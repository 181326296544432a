"""Per-cell semantics of computation strings on the GPU, in every kernel family: the programs of
``test_expr_lowering.py`` run on signed, seeded inputs with exact values planted at fixed cells.

Three tiers of reference:

* the table's compound strings against the oracle (``reference_numpy``), at the suite's tolerances;
* operations IEEE arithmetic rounds correctly (unary minus, fabs, min, max, floor, ceil, sqrt, the four
  arithmetic operators, selection, comparisons stored as 1.0 / 0.0): bit for bit against numpy in the field
  type, subnormal operands and results included -- a flush-to-zero or fast-math build fails here;
* transcendental functions: in ulps of the result, against numpy evaluated in float64 (float32 kernels) or in
  the 80-bit ``np.longdouble`` (float64 kernels) and rounded to the field type.

The cluster kernels share the one-operator kernels' cell code and must match them bit for bit."""
import json
import os
import zlib

import numpy as np
import pytest

import test_expr_lowering as tl

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-12}
# largest error in ulps each function may have: one above the maximum measured on a B200 (1000 W power limit;
# CUDA 12.9 NVRTC without fast math) over these inputs in every configuration, which was
# float32: sin 1, cos 1, tan 3, sinh 3, cosh 2, tanh 2, exp 2, log 1, pow 1, pow of negative bases 1;
# float64: sin 1, cos 1, tan 2, sinh 1, cosh 1, tanh 1, exp 1, log 1, pow 1, pow of negative bases 1
ULP_BOUND = {
    "float32": {"sin": 2, "cos": 2, "tan": 4, "sinh": 4, "cosh": 3, "tanh": 3, "exp": 3, "log": 2, "pow": 2,
                "powi": 2},
    "float64": {"sin": 2, "cos": 2, "tan": 3, "sinh": 2, "cosh": 2, "tanh": 2, "exp": 2, "log": 2, "pow": 2,
                "powi": 2},
}
TABLE_PROGRAMS = [n for n, (g, _) in tl.PROGRAMS.items() if g in tl.SCALAR]


@pytest.fixture(scope="module")
def gpu(native_lib):
    from stencilflow_b200 import runtime
    return runtime.Runtime.get()


def _planted(dt):
    """Integers, half-integers and their negatives, signed zeros, subnormals and the smallest normal."""
    fi = np.finfo(dt)
    sub, tiny = fi.smallest_subnormal, fi.tiny
    return np.array([0.0, -0.0, 0.5, -0.5, 1.0, -1.0, 1.5, -1.5, 2.0, -2.0, 0.25, -1.75, sub, -sub, 3 * sub, -3 * sub,
                     tiny / 2, -tiny / 4, tiny, -1.5 * tiny], dtype=dt)


def _plant(a, b, dt):
    """At runs of cells at the start, in the middle and at the end of the grid: ``a`` takes each planted value in
    two k-neighbouring cells; ``b`` equals ``a`` at the first (-a at the second, so sums and differences of
    subnormals are subnormal), except where that would divide zero by zero."""
    vals = _planted(dt)
    fa, fb = a.reshape(-1), b.reshape(-1)
    n = fa.size
    for base in (0, n // 3, 2 * n // 3, n - 3 * len(vals)):
        for q, v in enumerate(vals):
            c = base + 3 * q
            fa[c] = fa[c + 1] = v
            if fb is not None:
                fb[c], fb[c + 1] = (v, -v) if v != 0 else (dt(0.5), dt(-0.5))


def _positive(rng, shape, dt):
    p = rng.uniform(0.1, 4.0, size=shape).astype(dt)
    fi = np.finfo(dt)
    flat = p.reshape(-1)
    for q, v in enumerate((fi.smallest_subnormal, 3 * fi.smallest_subnormal, fi.tiny / 2, fi.tiny, 1.0, 4.0, 0.25)):
        flat[7 * q] = flat[flat.size // 2 + q] = v
    return p


def make_inputs(name, case):
    _, dtype, shape = case
    dt = np.dtype(dtype).type
    group = tl.PROGRAMS[name][0]
    # seeded by program, type and grid, not by configuration: the cluster run gets the one-operator run's inputs
    rng = np.random.default_rng(zlib.crc32("{}/{}/{}".format(name, dtype, shape).encode()))
    out = {}
    if group in ("signed", "exact"):
        out["a"] = rng.uniform(-2.0, 2.0, size=shape).astype(dt)
        out["b"] = rng.uniform(-2.0, 2.0, size=shape).astype(dt)
        _plant(out["a"], out["b"], dt)
    elif group == "positive":
        out["a"] = _positive(rng, shape, dt)
        out["b"] = _positive(rng, shape, dt)
    elif group == "pow":
        out["a"] = rng.uniform(0.5, 2.0, size=shape).astype(dt)              # bases (also of t)
        out["b"] = rng.integers(-3, 4, size=shape).astype(dt)                # integer exponents of negative bases
    if group == "exact":
        out["p"] = _positive(rng, shape, dt)
    if group == "transcendental":
        out["a"] = rng.uniform(-2.0, 2.0, size=shape).astype(dt)
        _plant(out["a"], np.zeros_like(out["a"]), dt)
        out["p"] = _positive(rng, shape, dt)
        out["q"] = rng.uniform(0.5, 2.0, size=shape).astype(dt)
        out["e"] = rng.uniform(-2.0, 2.0, size=shape).astype(dt)
        out["n"] = -rng.uniform(0.5, 2.0, size=shape).astype(dt)
        out["m"] = rng.integers(-3, 4, size=shape).astype(dt)
    if group in tl.SCALAR:
        out["s"] = dt(tl.SCALAR[group])
    return out


def _run(path, inputs, case, specialize=None):
    from oracle import reference_numpy as rn
    from stencilflow_b200.cuda_program import CudaProgram
    prog = CudaProgram(path, plan_options=tl.plan_options(case, path), specialize_scalars=specialize)
    try:
        tl.check_families(prog.plan, case)
        info = rn.ProgramInfo(rn.load_program(path))
        outs = {o: np.zeros(info.shape, dtype=info.field_type(o)) for o in info.outputs}
        args = {(k + "_host" if np.ndim(v) > 0 else k): v for k, v in inputs.items()}
        args.update({k + "_host": v for k, v in outs.items()})
        prog(**args)
    finally:
        prog.close()
    return outs


def _reference(path, inputs):
    from oracle import reference_numpy as rn
    with np.errstate(all="ignore"):
        return rn.run_reference(path, inputs)


def _trim(arr, halo):
    from oracle import reference_numpy as rn
    return rn.trim_halo(arr, halo)


def _run_case(name, case, tmp_path, monkeypatch, specialize=None):
    tl.clean_environment(monkeypatch, case)
    path, halos = tl.write_program(name, case, tmp_path)
    inputs = make_inputs(name, case)
    return path, halos, inputs, _run(path, inputs, case, specialize)


def _check_cluster_matches_general(name, case, tmp_path, monkeypatch, got, halos):
    if case[0] != "cluster":
        return
    general = ("general",) + tuple(case[1:])
    _, _, _, ref = _run_case(name, general, tmp_path, monkeypatch)
    for field, arr in got.items():
        assert _trim(arr, halos[field]).tobytes() == _trim(ref[field], halos[field]).tobytes(), field


def _check_oracle(path, halos, inputs, got, case):
    """At the suite's tolerances.  Inputs and results are of order one and cross zero, so near zero the bound is
    absolute at that scale: |got - ref| <= tol * max(|ref|, 1)."""
    expected = _reference(path, inputs)
    for field, ref in expected.items():
        r = _trim(ref, halos[field]).astype(np.float64)
        g = _trim(got[field], halos[field]).astype(np.float64)
        assert np.isfinite(r).all(), field
        err = np.abs(r - g) / np.maximum(np.abs(r), 1.0)
        worst = np.unravel_index(np.nanargmax(np.where(np.isnan(err), np.inf, err)), err.shape)
        assert np.isfinite(g).all() and err.max() <= TOL[case[1]], \
            "{} {}: err {} at {}: got {} want {}".format(tl.case_id(case), field, err[worst], worst, g[worst], r[worst])


@pytest.mark.parametrize("name", TABLE_PROGRAMS)
@pytest.mark.parametrize("case", tl.CASES, ids=tl.case_id)
def test_table_matches_the_oracle(gpu, tmp_path, monkeypatch, case, name):
    path, halos, inputs, got = _run_case(name, case, tmp_path, monkeypatch)
    _check_oracle(path, halos, inputs, got, case)
    _check_cluster_matches_general(name, case, tmp_path, monkeypatch, got, halos)


@pytest.mark.parametrize("name", TABLE_PROGRAMS)
@pytest.mark.parametrize("case", [c for c in tl.CASES if c[2] == tl.SMALL and c[0] in ("general", "packed", "stream64")],
                         ids=tl.case_id)
def test_specialized_scalars_match_the_oracle(gpu, tmp_path, monkeypatch, case, name):
    """``s`` as a literal of the kernel (the compiler may then fold and contract differently, so not bit for bit
    the kernel with ``s`` as a parameter)."""
    group = tl.PROGRAMS[name][0]
    path, halos, inputs, got = _run_case(name, case, tmp_path, monkeypatch, specialize={"s": tl.SCALAR[group]})
    _check_oracle(path, halos, inputs, got, case)


@pytest.mark.parametrize("case", tl.CASES, ids=tl.case_id)
def test_correctly_rounded_operations_are_exact(gpu, tmp_path, monkeypatch, case):
    path, halos, inputs, got = _run_case("exact", case, tmp_path, monkeypatch)
    dt = np.dtype(case[1]).type
    # numpy in the field type, with subnormals (copy boundaries keep the oracle there)
    expected = _reference(path, inputs)
    fi = np.finfo(dt)
    a = inputs["a"]
    assert ((np.abs(a) < fi.tiny) & (a != 0)).sum() >= 16
    bad = []
    for field, ref in expected.items():
        assert ref.dtype == dt
        if not np.array_equal(ref, got[field]):
            diff = np.argwhere(ref != got[field])
            c = tuple(diff[0])
            bad.append("{}: {} cells, first {} got {!r} want {!r}".format(field, len(diff), c, got[field][c], ref[c]))
    # subnormal results survive
    sub = (np.abs(expected["min"]) < fi.tiny) & (expected["min"] != 0)
    assert sub.any()
    assert not bad, bad
    _check_cluster_matches_general("exact", case, tmp_path, monkeypatch, got, halos)


def _ulps(got, ref):
    """|got - ref| in units of the last place of ``ref`` (both of the field type)."""
    ref64 = ref.astype(np.float64)
    return np.abs(got.astype(np.float64) - ref64) / np.spacing(np.abs(ref)).astype(np.float64)


def test_ulps_of_correctly_rounded_values():
    x = np.float32(1.5)
    assert _ulps(np.array([np.nextafter(x, np.float32(2))]), np.array([x]))[0] == 1.0
    sub = np.finfo(np.float64).smallest_subnormal
    assert _ulps(np.array([3 * sub]), np.array([sub]))[0] == 2.0


@pytest.mark.parametrize("case", tl.CASES, ids=tl.case_id)
def test_transcendental_functions_within_their_ulp_bounds(gpu, tmp_path, monkeypatch, case):
    path, halos, inputs, got = _run_case("transcendental", case, tmp_path, monkeypatch)
    dtype = case[1]
    dt = np.dtype(dtype).type
    wide = np.float64 if dtype == "float32" else np.longdouble
    x = {k: v.astype(wide) for k, v in inputs.items()}
    exact = {"sin": np.sin(x["a"]), "cos": np.cos(x["a"]), "tan": np.tan(x["a"]), "sinh": np.sinh(x["a"]),
             "cosh": np.cosh(x["a"]), "tanh": np.tanh(x["a"]), "exp": np.exp(x["a"]), "log": np.log(x["p"]),
             "pow": np.power(x["q"], x["e"]), "powi": np.power(x["n"], x["m"])}
    measured, bad = {}, []
    for fn, want in exact.items():
        ref = want.astype(dt)
        assert np.isfinite(ref).all() and np.isfinite(got[fn]).all(), fn
        ulps = _ulps(got[fn], ref)
        measured[fn] = float(ulps.max())
        if measured[fn] > ULP_BOUND[dtype][fn]:
            c = np.unravel_index(np.argmax(ulps), ulps.shape)
            bad.append("{}: {} ulp at {}: x={!r} got {!r} want {!r}".format(fn, measured[fn], c,
                                                                         [inputs[k][c] for k in ("a", "p", "q", "e", "n", "m")],
                                                                         got[fn][c], ref[c]))
    print("ulp maxima", tl.case_id(case), measured)
    assert not bad, bad
    _check_cluster_matches_general("transcendental", case, tmp_path, monkeypatch, got, halos)


@pytest.mark.parametrize("unroll", ["1", "6"])
def test_copy_boundaries_on_a_grid_with_boundary_free_trips(gpu, tmp_path, monkeypatch, unroll):
    """The copy-boundary Jacobi-3D chain of the test programs on a grid whose fused pass runs trips without boundary
    code: the last operator's i-1 tap at plane 0 must read its own plane, not one outside the domain.  Against the
    oracle and, bit for bit, the one-operator kernels."""
    from conftest import program_path
    from oracle import reference_numpy as rn
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    for k in [k for k in os.environ if k.startswith("SFB200_") and k != "SFB200_CACHE"]:
        monkeypatch.delenv(k)
    monkeypatch.setenv("SFB200_UNROLL", unroll)
    with open(program_path("jacobi3d_12x12x16_3itr_copy")) as f:
        desc = json.load(f)
    shape = [24, 200, 384]
    desc["dimensions"] = shape
    path = str(tmp_path / "jacobi3d_copy_large.json")
    with open(path, "w") as f:
        json.dump(desc, f)
    a = np.random.default_rng(3).uniform(0.0, 1.0, size=shape).astype(np.float32)
    expected = rn.run_reference(path, {"a": a})["b2"]
    results = {}
    for label, opts in (("unfused", PlanOptions(fuse=False)), ("fused", PlanOptions(max_depth=3))):
        prog = CudaProgram(path, plan_options=opts)
        try:
            streamed = [l for l in prog.lowered.launches if l.family == "streamed"]
            if label == "fused":
                assert len(streamed) == 1
                rows, cols = streamed[0].info["tile"]
                assert shape[1] >= 3 * rows and shape[2] >= 3 * cols
            out = np.zeros(shape, np.float32)
            prog(a_host=a, b2_host=out)
        finally:
            prog.close()
        err = rn.max_relative_error(expected, out)
        assert err <= TOL["float32"], "{}: max rel err {} at {}".format(
            label, err, np.unravel_index(np.argmax(np.abs(expected - out)), shape))
        results[label] = out.tobytes()
    assert results["fused"] == results["unfused"]

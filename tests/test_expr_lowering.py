"""Computation strings through every per-cell emitter (no GPU): a table of strings that covers the grammar of
``expr.py``, lowered in each kernel family and compiled with NVRTC.  ``test_expr_semantics_gpu.py`` runs the same
programs on the GPU against the oracle.

Each table string is the consumer of an intermediate ``t = a[i,j,k]``, so that in a fused pass it reads ``t``
through the exchange ring; its taps reach the i, j and k boundaries under constant, shrink and copy conditions.
Independent consumers of one producer share a program to keep the number of compiles down."""
import json
import os
import re

import pytest


DIMS = ["i", "j", "k"]
SCALAR = {"signed": -0.75, "positive": 1.25, "pow": 1.5}     # the 0-D input ``s`` of each input group
C0 = 0.25                                                     # the program constant ``c0``

# (consumer name, input group, computation string).  The groups fix the input ranges (test_expr_semantics_gpu):
# "signed" [-2, 2], "positive" [0.1, 4] (log, sqrt), "pow" bases in [0.5, 2] and integer-valued exponents.
# Literals the float32 and float64 lowerings could round differently are kept dyadic.
TABLE = [
    ("trig", "signed",
     "r = sin(t[i-1,j,k]) + cos(t[i,j+1,k]) * tan(0.5 * a[i,j,k-1]) - sin(s) * cos(t[i,j,k])"),
    ("hyper", "signed",
     "r = sinh(t[i,j,k]) - cosh(a[i+1,j,k]) * 0.25 + tanh(t[i,j-1,k+1] * s) + tanh(c0)"),
    ("expround", "signed",
     "r = exp(t[i,j,k-1]) * 0.25 + floor(t[i+1,j,k] * 4.0) - ceil(b[i,j+1,k] * 2.0) + floor(t[i,j,k]) "
     "+ ceil(a[i,j,k]) + fabs(t[i,j,k+1]) - abs(a[i,j,k]) + abs(s) + exp(c0)"),
    ("minmax", "signed",
     "r = min(t[i,j,k], s) + max(c0, a[i,j+1,k]) + min(a[i-1,j,k], t[i,j,k+1]) + max(t[i,j,k-1], b[i,j,k]) "
     "+ min(s, c0) + max(b[i,j,k], s)"),
    ("compare", "signed",
     "r = (1.0 if t[i,j,k] < a[i,j,k+1] else 0.0) + (2.0 if t[i-1,j,k] <= 0.5 else 0.0) "
     "+ (4.0 if t[i,j+1,k] > b[i,j,k] else 0.0) + (8.0 if a[i,j,k+1] >= -0.25 else 0.0) "
     "+ (16.0 if t[i,j,k] == b[i,j,k] else 0.0) + (32.0 if t[i,j,k-1] != a[i,j,k] else 0.0) "
     "+ (64.0 if s < c0 else 0.0)"),
    ("logic", "signed",
     "c = t[i,j,k] > 0.5 and a[i,j-1,k] < 0.25 and b[i,j,k] > -0.5; "
     "d = t[i+1,j,k] < -0.5 or a[i,j,k] > 1.5 or not (b[i,j,k+1] <= 0.25); "
     "e = not (s > c0) or t[i,j,k] == a[i,j,k]; "
     "r = (1.0 if c else 0.0) + (2.0 if d else 0.0) + (4.0 if not c else 0.0) + (8.0 if e else 0.0)"),
    ("select", "signed",
     "c = (t[i,j,k] > 0.5) if a[i,j,k] > 0.0 else (t[i,j,k-1] < 0.25); "
     "r = t[i,j,k] if c else (b[i-1,j,k] if t[i,j+1,k] < 0.0 else (-a[i,j,k] if s > c0 else 2.0))"),
    ("negate", "signed",
     "x = t[i,j,k] * 0.5; y = -s; r = -t[i-1,j,k] + y * a[i,j,k-1] - (-x) + -(c0 * s) - -b[i,j+1,k]"),
    # the FMA shapes of the packed emitter, the uniform operand in each position it can take; the odd k-offsets
    # are not register pairs and take the conventional path
    ("fma_add", "signed",
     "p1 = s * t[i,j,k] + a[i,j,k]; p2 = t[i,j,k] * s + b[i,j,k]; p3 = t[i,j,k] * a[i,j,k] + c0; "
     "p4 = t[i,j,k] * a[i,j,k] + b[i,j,k]; p5 = a[i,j,k] + s * t[i,j,k]; p6 = b[i,j,k] + t[i,j,k] * c0; "
     "p7 = s + t[i,j,k] * b[i,j,k]; p8 = t[i-1,j,k] + t[i,j,k+1] * a[i,j+1,k]; "
     "r = p1 + p2 + p3 + p4 + p5 + p6 + p7 + p8"),
    ("fma_sub", "signed",
     "m1 = t[i,j,k] * a[i,j,k] - s; m2 = s * t[i,j,k] - b[i,j,k]; m3 = t[i,j,k] * c0 - a[i,j,k]; "
     "m4 = t[i,j,k] * a[i,j,k] - b[i,j-1,k]; n1 = s - t[i,j,k] * b[i,j,k]; n2 = a[i,j,k] - c0 * t[i,j,k]; "
     "n3 = b[i,j,k] - t[i,j,k] * s; n4 = b[i+1,j,k] - t[i,j,k] * a[i,j,k-1]; "
     "r = m1 + 2.0 * m2 + 4.0 * m3 + 8.0 * m4 + 0.5 * n1 + 0.25 * n2 - n3 - 2.0 * n4"),
    ("uniform_temps", "signed",
     "u = s * c0; v = u + 2.0; w = -u; z = 3.0; "
     "r = t[i,j,k] * v + (u if s > c0 else w) + a[i,j+1,k] * w - z * t[i,j,k-1] + b[i-1,j,k]"),
    ("reassign", "signed",
     "x = t[i,j,k]; x = x + t[i,j,k+1]; x = x * 0.5; y = a[i-1,j,k]; y = y - x; r = x - y * b[i,j+1,k]"),
    ("bool_reassign", "signed",
     "c = t[i,j,k] > 0.5; c = c and a[i,j,k] < 0.75; c = c or b[i,j+1,k] < -1.5; "
     "r = 1.0 if c else 2.0 + t[i-1,j,k-1]"),
    ("retype", "signed",
     "c = t[i,j,k] > 0.5; c = t[i,j,k] * 2.0 + a[i+1,j,k]; d = t[i,j,k] * 2.0; d = d > a[i,j-1,k]; "
     "r = c + d + (1.0 if d else -1.0) - t[i,j,k+1]"),
    # the result is the last statement's target, not the operator's name
    ("named", "signed",
     "x = t[i,j,k] + a[i,j,k+1]; y = x * x - b[i-1,j,k] + t[i,j-1,k]"),
    ("literals", "signed",
     "r = t[i,j,k] * 1e-3 + 2 * a[i,j,k] + (1 / 2) * b[i,j-1,k] + (1.0 if True else 0.0) + 3 "
     "+ (0.5 if False else t[i+1,j,k]) - 1.5e1 * c0 + t[i,j,k+1]"),
    ("logsqrt", "positive",
     "r = log(t[i,j,k]) + sqrt(a[i,j+1,k]) * log(b[i-1,j,k]) - sqrt(t[i,j,k-1] * s) + log(s) + sqrt(c0)"),
    ("powers", "pow",
     "r = pow(t[i,j,k], s) + pow(a[i,j+1,k], t[i,j,k-1]) + pow(-t[i-1,j,k], 3.0) + pow(-t[i,j,k], b[i,j,k]) "
     "+ pow(c0, t[i,j,k+1]) + pow(s, c0)"),
]

# operations that are correctly rounded in IEEE arithmetic: one operator each, no literal, copy boundaries only
# (they keep the oracle in the field type), compared bit for bit
EXACT = [
    ("neg", "-a[i,j,k]"), ("fabs", "fabs(a[i,j,k])"), ("abs", "abs(b[i,j,k])"),
    ("min", "min(a[i,j,k], b[i,j,k])"), ("max", "max(a[i,j,k], b[i,j,k])"),
    ("floor", "floor(a[i,j,k])"), ("ceil", "ceil(b[i,j,k])"), ("sqrt", "sqrt(p[i,j,k])"),
    ("add", "a[i,j,k] + b[i,j,k]"), ("sub", "a[i,j,k] - b[i,j,k]"), ("mul", "a[i,j,k] * b[i,j,k]"),
    ("div", "a[i,j,k] / b[i,j,k]"), ("subk", "a[i,j,k+1] - a[i,j,k]"), ("addj", "b[i,j-1,k] + b[i,j,k]"),
    ("sel", "a[i,j,k] if a[i,j,k] < b[i,j,k] else b[i,j,k]"),
    ("lt", "a[i,j,k] < b[i,j,k]"), ("le", "a[i,j,k] <= b[i,j,k]"), ("gt", "a[i,j,k] > b[i,j,k]"),
    ("ge", "a[i,j,k] >= b[i,j,k]"), ("eq", "a[i,j,k] == b[i,j,k]"), ("ne", "a[i,j,k] != b[i,j,k]"),
]

# transcendental functions, one operator each, measured in ulps of the result
TRANSCENDENTAL = [
    ("sin", "sin(a[i,j,k])"), ("cos", "cos(a[i,j,k])"), ("tan", "tan(a[i,j,k])"), ("sinh", "sinh(a[i,j,k])"),
    ("cosh", "cosh(a[i,j,k])"), ("tanh", "tanh(a[i,j,k])"), ("exp", "exp(a[i,j,k])"), ("log", "log(p[i,j,k])"),
    ("pow", "pow(q[i,j,k], e[i,j,k])"), ("powi", "pow(n[i,j,k], m[i,j,k])"),
]

SMALL = [12, 20, 32]
# float32 / float64 grids on which the fused passes have tiles whose halo lies inside the domain (boundary-free trips)
LARGE = {"float32": [20, 200, 384], "float64": [20, 200, 256]}
UNALIGNED = {"float32": [12, 20, 30], "float64": [12, 20, 31]}   # innermost rows of 120 and 248 bytes

# label -> (PlanOptions keywords, environment, intended family); max_depth None = as many as the program has.
# The fused passes are not unrolled over streamed steps: the cell code is the same, the source a sixth as long
# (NVRTC time dominates these tests).
ONE_STEP = {"SFB200_UNROLL": "1"}
CONFIGS = {
    "general": (dict(fuse=False), {}, "general"),
    "packed": (dict(max_depth=None), ONE_STEP, "streamed"),
    "scalar": (dict(max_depth=None), dict(ONE_STEP, SFB200_PACK="0"), "streamed"),
    "stream64": (dict(max_depth=None), ONE_STEP, "streamed"),
    "unaligned": (dict(max_depth=None, unaligned=1), ONE_STEP, "streamed"),
    "cluster": (dict(cluster=1), {}, "cluster"),
}
# (configuration, dtype, shape)
CASES = [
    ("general", "float32", SMALL), ("general", "float64", SMALL),
    ("packed", "float32", SMALL), ("packed", "float32", LARGE["float32"]),
    ("scalar", "float32", SMALL),
    ("stream64", "float64", SMALL), ("stream64", "float64", LARGE["float64"]),
    ("unaligned", "float32", UNALIGNED["float32"]), ("unaligned", "float64", UNALIGNED["float64"]),
    ("cluster", "float32", SMALL), ("cluster", "float64", SMALL),
]
CONSUMERS_PER_PROGRAM = 5


def case_id(case):
    config, dtype, shape = case
    return "{}-{}-{}".format(config, dtype, "x".join(map(str, shape)))


def _groups():
    """Table programs: (name, group, [(consumer, string)]), at most CONSUMERS_PER_PROGRAM consumers each."""
    out = []
    for group in SCALAR:
        rows = [(n, cs) for n, g, cs in TABLE if g == group]
        for p in range(0, len(rows), CONSUMERS_PER_PROGRAM):
            out.append(("{}{}".format(group, p // CONSUMERS_PER_PROGRAM), group, rows[p:p + CONSUMERS_PER_PROGRAM]))
    return out


PROGRAMS = {name: (group, rows) for name, group, rows in _groups()}
PROGRAMS["exact"] = ("exact", [(n, "{} = {}".format(n, cs)) for n, cs in EXACT])
PROGRAMS["transcendental"] = ("transcendental", [(n, "{} = {}".format(n, cs)) for n, cs in TRANSCENDENTAL])

INPUTS = {"signed": ["a", "b"], "positive": ["a", "b"], "pow": ["a", "b"],
          "exact": ["a", "b", "p"], "transcendental": ["a", "p", "q", "e", "n", "m"]}


def parse(cs):
    from stencilflow_b200 import expr
    dims = {f: list(DIMS) for f in ("t", "a", "b", "p", "q", "e", "n", "m")}
    dims["s"] = []
    return expr.parse_computation(cs, dims, DIMS)


def _boundaries(cs, n):
    """Boundary conditions of consumer ``n``: constant, shrink and copy rotate over t, a and b (copy only where
    the centre tap is read, which a copy boundary needs).  Returns (conditions, halo to trim)."""
    from stencilflow_b200 import expr
    kinds = ("constant", "shrink", "copy")
    taps = expr.collect_taps(parse(cs))
    bcs, halo = {}, 0
    for m, field in enumerate(sorted(taps)):
        offsets = taps[field]
        if not any(any(o) for o in offsets):
            continue
        kind = kinds[(n + m) % 3]
        if kind == "copy" and (0, 0, 0) not in offsets:
            kind = "constant"
        bcs[field] = {"type": "copy"} if kind == "copy" else (
            {"type": "shrink"} if kind == "shrink" else {"type": "constant", "value": 0.5})
        if kind == "shrink":
            halo = max([halo] + [abs(o) for off in offsets for o in off])
    return bcs, halo


def program_desc(name, dtype, shape):
    """JSON description of table program ``name`` and {output: halo}."""
    from stencilflow_b200 import expr
    group, rows = PROGRAMS[name]
    inputs = {f: {"data": "constant:0.5", "data_type": dtype} for f in INPUTS[group]}
    ops, halos = {}, {}
    if group in SCALAR:
        inputs["s"] = {"data": SCALAR[group], "data_type": dtype, "input_dims": []}
        ops["t"] = {"computation_string": "t = a[i,j,k]", "data_type": dtype, "boundary_conditions": {}}
        for n, (consumer, cs) in enumerate(rows):
            bcs, halos[consumer] = _boundaries(cs, n)
            ops[consumer] = {"computation_string": cs, "data_type": dtype, "boundary_conditions": bcs}
    else:
        for consumer, cs in rows:
            fields = {f for f, offs in expr.collect_taps(parse(cs)).items() if any(any(o) for o in offs)}
            ops[consumer] = {"computation_string": cs, "data_type": dtype,
                             "boundary_conditions": {f: {"type": "copy"} for f in sorted(fields)}}
            halos[consumer] = 0
    desc = {"inputs": inputs, "outputs": [o for o in ops if o != "t"], "dimensions": list(shape), "program": ops}
    if group in SCALAR:
        desc["constants"] = {"c0": {"data_type": dtype, "value": C0}}
    return desc, halos


def write_program(name, case, directory):
    config, dtype, shape = case
    desc, halos = program_desc(name, dtype, shape)
    path = os.path.join(str(directory), "{}_{}.json".format(name, case_id(case)))
    with open(path, "w") as f:
        json.dump(desc, f)
    return path, halos


def plan_options(case, path):
    from stencilflow_b200.planner import PlanOptions
    opts = dict(CONFIGS[case[0]][0])
    if "max_depth" in opts:
        with open(path) as f:
            opts["max_depth"] = len(json.load(f)["program"])
    return PlanOptions(**opts)


def clean_environment(monkeypatch, case):
    for k in list(os.environ):
        if k.startswith("SFB200_") and k != "SFB200_CACHE":
            monkeypatch.delenv(k)
    for k, v in CONFIGS[case[0]][1].items():
        monkeypatch.setenv(k, v)


def check_families(plan, case):
    """The launches are of the family the configuration is for."""
    config, dtype, shape = case
    family = CONFIGS[config][2]
    launches = plan.lowered.launches
    assert launches and all(l.family == family for l in launches), [l.family for l in launches]
    if family == "cluster":
        assert len(launches) == 1
    if config == "unaligned":
        assert all(l.info.get("unaligned") for l in launches)
    if shape == LARGE.get(dtype) and family == "streamed":
        for l in launches:
            rows, cols = l.info["tile"]
            assert shape[1] >= 3 * rows and shape[2] >= 3 * cols, (l.info["tile"], shape)


def _lower(name, case, tmp_path, monkeypatch, specialize=None):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.planner import plan_program
    from stencilflow_b200.stencil_op import make_program
    clean_environment(monkeypatch, case)
    path, _ = write_program(name, case, tmp_path)
    plan = plan_program(make_program(KernelChainGraph(path)), plan_options(case, path), specialize=specialize)
    check_families(plan, case)
    return path, plan


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_table_lowers_to_the_family_and_compiles(native_lib, tmp_path, monkeypatch, case):
    from stencilflow_b200.cuda_program import CudaProgram
    monkeypatch.setenv("SFB200_CACHE", str(tmp_path / "cache"))
    for name in PROGRAMS:
        path, plan = _lower(name, case, tmp_path, monkeypatch)
        prog = CudaProgram(path, plan_options=plan_options(case, path), allocate=False)
        assert len(prog.image) > 0, name
        assert prog.lowered.source == plan.lowered.source, name


@pytest.mark.parametrize("case", [c for c in CASES if c[2] == SMALL and c[0] in ("general", "packed", "stream64")],
                         ids=case_id)
def test_specialized_scalars_compile(native_lib, tmp_path, monkeypatch, case):
    """The 0-D input as a literal of the kernel (``specialize_scalars``) rather than a kernel parameter."""
    from stencilflow_b200.cuda_program import CudaProgram
    monkeypatch.setenv("SFB200_CACHE", str(tmp_path / "cache"))
    for name, (group, _) in PROGRAMS.items():
        if group not in SCALAR:
            continue
        path, plan = _lower(name, case, tmp_path, monkeypatch, specialize={"s": SCALAR[group]})
        assert not [a for l in plan.lowered.launches for a in l.args if a[0] == "scalar"], name
        prog = CudaProgram(path, plan_options=plan_options(case, path), specialize_scalars={"s": SCALAR[group]},
                           allocate=False)
        assert len(prog.image) > 0, name


@pytest.mark.parametrize("string", [
    "c = t[i,j,k] > 0.5; c = c and a[i,j,k] < 0.7; r = 1.0 if c else 2.0",
    "x = t[i,j,k]; x = x + t[i,j,k+1]; x = x * 0.5; r = x",
])
@pytest.mark.parametrize("case", [c for c in CASES if c[2] == SMALL or c[0] == "unaligned"], ids=case_id)
def test_reassigned_temporaries_compile(native_lib, tmp_path, monkeypatch, case, string):
    """Two strings that once failed to compile: a boolean temporary assigned twice (an assignment to a const
    bool) in the one-operator and cluster kernels, and a temporary assigned three times (a name declared
    twice) in the float64 and one-cell-at-a-time fused passes."""
    from stencilflow_b200.cuda_program import CudaProgram
    monkeypatch.setenv("SFB200_CACHE", str(tmp_path / "cache"))
    clean_environment(monkeypatch, case)
    config, dtype, shape = case
    desc = {"inputs": {"a": {"data": "constant:0.5", "data_type": dtype}}, "outputs": ["r"],
            "dimensions": list(shape),
            "program": {"t": {"computation_string": "t = a[i,j,k]", "data_type": dtype, "boundary_conditions": {}},
                        "r": {"computation_string": string, "data_type": dtype,
                              "boundary_conditions": {"t": {"type": "constant", "value": 0.0}}}}}
    path = str(tmp_path / "reassign.json")
    with open(path, "w") as f:
        json.dump(desc, f)
    prog = CudaProgram(path, plan_options=plan_options(case, path), allocate=False)
    check_families(prog.plan, case)
    assert len(prog.image) > 0


def test_reassignment_takes_the_type_of_its_own_value():
    """A number assigned to a name that held a boolean stays a number (and the reverse), in every emitter that
    declares C variables."""
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.planner import PlanOptions, plan_program
    from stencilflow_b200.stencil_op import make_program
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        path, _ = write_program("signed2", ("general", "float64", SMALL), d)
        src = plan_program(make_program(KernelChainGraph(path)), PlanOptions(fuse=False)).lowered.source
    # retype: c bool then double, d double then bool
    assert re.search(r"const bool v0_t(\d+) = .*\n  double v0_t\1_1 = ", src)
    assert re.search(r"  double v0_t(\d+) = .*\n(  .*\n)*?  const bool v0_t\1_1 = ", src)


def _constructs(stmts):
    from stencilflow_b200 import expr as ex
    seen = set()
    for s in stmts:
        for e in ex.walk(s.value):
            if isinstance(e, ex.Call):
                seen.add(("call", e.fn))
                if len(e.args) == 2:
                    kinds = {"field" if any(isinstance(x, ex.Tap) for x in ex.walk(a)) else "uniform" for a in e.args}
                    if kinds == {"field", "uniform"}:
                        seen.add(("mixed call", e.fn))
            elif isinstance(e, ex.Cmp):
                seen.add(("cmp", e.op))
            elif isinstance(e, ex.Logic):
                seen.add(("logic", e.op, min(len(e.args), 3)))
            elif isinstance(e, ex.Select):
                seen.add("select")
                if isinstance(e.a, ex.Select) or isinstance(e.b, ex.Select):
                    seen.add("nested select")
                if all(isinstance(x, (ex.Cmp, ex.Logic)) for x in (e.a, e.b)):
                    seen.add("boolean select")
            elif isinstance(e, ex.Neg):
                seen.add(("neg", type(e.a).__name__))
            elif isinstance(e, ex.Const):
                seen.add(("literal", type(e.value).__name__))
    return seen


def test_table_covers_the_grammar():
    """Every function (both spellings of fabs), comparison, logic operator, ternary shape and literal kind appears
    in the table: a function or operator added to ``expr.py`` without a case here fails this test."""
    from stencilflow_b200 import expr as ex
    seen = set()
    for _, _, cs in TABLE:
        seen |= _constructs(parse(cs))
    need = {("call", f) for f in ex.FUNCTIONS}
    need |= {("mixed call", f) for f, (_, arity) in ex.FUNCTIONS.items() if arity == 2}
    need |= {("cmp", op) for op in ex._CMPOPS.values()}
    need |= {("logic", "and", 3), ("logic", "or", 3), ("logic", "not", 1)}
    need |= {"select", "nested select", "boolean select"}
    need |= {("neg", "Tap"), ("neg", "Var"), ("neg", "Bin")}
    need |= {("literal", "int"), ("literal", "float"), ("literal", "bool")}
    assert need <= seen, sorted(map(str, need - seen))
    strings = [cs for _, _, cs in TABLE]
    assert any("1e-3" in cs for cs in strings) and any("(1 / 2)" in cs for cs in strings)
    # the exact and transcendental programs cover their functions too
    exact = set().union(*(_constructs(parse("r = " + cs)) for _, cs in EXACT))
    assert {("call", f) for f in ("fabs", "abs", "min", "max", "floor", "ceil", "sqrt")} <= exact
    assert {("cmp", op) for op in ex._CMPOPS.values()} <= exact
    trans = set().union(*(_constructs(parse("r = " + cs)) for _, cs in TRANSCENDENTAL))
    assert {("call", f) for f in ("sin", "cos", "tan", "sinh", "cosh", "tanh", "exp", "log", "pow")} <= trans


def test_table_temporaries():
    """Temporaries from uniform values only, assigned two and three times, booleans reassigned, reassignments that
    change the type both ways, and a result named other than its operator."""
    stmts = {n: parse(cs) for n, _, cs in TABLE}
    counts = {n: {t: [s.target for s in st].count(t) for t in {s.target for s in st}} for n, st in stmts.items()}
    assert any(3 in c.values() for c in counts.values()) and any(2 in c.values() for c in counts.values())
    from stencilflow_b200 import expr as ex

    def is_bool(e):
        return isinstance(e, (ex.Cmp, ex.Logic))
    changes = set()
    for st in stmts.values():
        last = {}
        for s in st:
            if s.target in last:
                changes.add((last[s.target], is_bool(s.value)))
            last[s.target] = is_bool(s.value)
    assert {(True, True), (True, False), (False, True), (False, False)} <= changes
    assert any(not any(isinstance(e, ex.Tap) for e in ex.walk(s.value)) and
               any(isinstance(e, ex.Var) for e in ex.walk(s.value)) for st in stmts.values() for s in st)
    assert any(st[-1].target not in ("r",) for st in stmts.values())


def test_every_consumer_reaches_the_boundaries_under_each_condition():
    kinds = set()
    for name, (group, rows) in PROGRAMS.items():
        if group not in SCALAR:
            continue
        desc, _ = program_desc(name, "float32", SMALL)
        for consumer, cs in rows:
            from stencilflow_b200 import expr
            taps = expr.collect_taps(parse(cs))
            assert "t" in taps, consumer
            reach = [any(off[d] for offs in taps.values() for off in offs) for d in range(3)]
            assert all(reach), (consumer, reach)
            kinds |= {bc["type"] for bc in desc["program"][consumer]["boundary_conditions"].values()}
    assert kinds == {"constant", "shrink", "copy"}


def test_packed_emitter_branches(tmp_path, monkeypatch):
    """The float32 fused passes of the table together use every kind of value of the packed emitter: packed FMA,
    addition, subtraction and multiplication, a uniform operand widened to a pair, and boolean lane pairs."""
    sources = []
    for case in CASES:
        if case[0] != "packed":
            continue
        for name in PROGRAMS:
            sources.append(_lower(name, case, tmp_path, monkeypatch)[1].lowered.source)
    text = "\n".join(sources)
    for fn in ("sf_fma2(", "sf_add2(", "sf_sub2(", "sf_mul2("):
        assert fn in text, fn
    assert re.search(r"make_float2\(([^,]+), \1\)", text)
    assert re.search(r"const bool (\w+)l = \(.*\), \1h = \(", text)

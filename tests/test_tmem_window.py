"""Tensor-memory window slots of the fused 3-D pass (no GPU): which slots qualify, what the register estimate
and the shared-memory budget make of them, and what the generator emits."""
import pytest

from conftest import program_path


def _program(name):
    return _program_at(program_path(name))


def _program_at(path):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    return make_program(KernelChainGraph(path))


def _analysis(prog, ops=None):
    from stencilflow_b200 import lower_stream
    return lower_stream.GroupAnalysis(prog, ops or list(prog.ops), exchange_cols=False)


def _config1():
    from stencilflow_b200 import programs
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    name, prog, _ = programs.baseline_config(1)
    return make_program(KernelChainGraph(programs.write_program(prog, name)))


def test_jacobi3d_parks_the_oldest_plane_of_every_window():
    """A 7-point chain reads the i-1 plane of each window only at the consumer's own cell: all four windows
    of a 4-operator pass qualify, at age 2; the last result is not consumed and has no window."""
    prog = _program("ref_jacobi3d_32x32x32_8itr")
    ana = _analysis(prog, list(prog.ops)[:4])
    assert {n: i.window for n, i in ana.fields.items() if i.consumed} == {n: 3 for n in ana.tmem_ages}
    assert len(ana.tmem_ages) == 4 and set(ana.tmem_ages.values()) == {2}


def test_hdiff_parks_only_the_planes_read_at_the_own_cell():
    """hdiff streamed along i: the i+1 tap of ``lap`` makes ``inp`` four planes deep and ``flx`` three; their
    oldest planes are read at the own cell only.  ``lap`` and ``fly`` end on planes read by j-neighbours."""
    ana = _analysis(_program("hdiff_24x28x16"))
    assert dict(ana.tmem_ages) == {"inp": 3, "flx": 2}
    assert ana.fields["lap"].window == 2 and ana.fields["fly"].window == 2


@pytest.mark.parametrize("name", ["jacobi2d_64x64_4itr_const_f32", "jacobi2d_96x128_6itr_shrink_f64"])
def test_no_tensor_memory_in_2d_passes(name):
    """2-D passes run several CTAs per SM: whatever their windows, they never get tensor memory."""
    from stencilflow_b200 import lower_stream
    ana = _analysis(_program(name))
    built = 0
    for V in (2, 4):
        for (R, WR, WC, KS) in [(1, 1, 1, 32), (1, 1, 2, 32), (1, 1, 8, 32)]:
            try:
                geo = lower_stream.Geometry(ana, V, R, WR, WC, 2, KS, tmem=True)
            except lower_stream.NotStreamable:
                continue
            built += 1
            assert not geo.tmem and geo.tmem_cols == 0
    assert built


def test_register_estimate_drops_by_the_parked_planes():
    prog = _config1()
    ana = _analysis(prog, list(prog.ops)[:4])
    assert ana.register_estimate(3, 4) == 168
    assert ana.register_estimate(3, 4, tmem=True) == 168 - 4 * 12
    assert ana.register_estimate(4, 4, tmem=True) == ana.register_estimate(4, 4) - 4 * 16


def test_r4_geometry_fits_shared_memory_and_tensor_memory():
    """R = 4 x 12 warps (24 row groups of 16 threads, a 96 x 64 tile), TMA ring 4 ahead: 221 KB of shared memory,
    and registers only with the planes parked; 16-word planes, two per field, four fields = the 128 columns
    of each warp."""
    from stencilflow_b200 import lower_stream
    prog = _config1()
    ana = _analysis(prog, list(prog.ops)[:4])
    geo = lower_stream.Geometry(ana, 4, 4, 24, 1, 4, 16, tmem=True)
    assert geo.tmem and geo.tmem_cols == 16 and 2 * geo.tmem_cols * len(ana.tmem_ages) == 128
    assert geo.smem == 221320 <= lower_stream.SMEM_LIMIT
    assert lower_stream.resident_estimate(geo) == 1
    assert ana.register_estimate(4, 4, tmem=True) <= lower_stream.register_limit(geo.NT) < ana.register_estimate(4, 4)
    assert lower_stream.Geometry(ana, 4, 4, 24, 1, 4, 16).smem == geo.smem - 16


def test_generated_pass_allocates_parks_fetches_and_frees():
    from stencilflow_b200 import lower_stream
    prog = _config1()
    ops = list(prog.ops)[:4]
    ana = _analysis(prog, ops)
    geo = lower_stream.Geometry(ana, 4, 3, 24, 1, 5, 16, tmem=True)
    gen = lower_stream.StreamKernelGen(prog, ops, ana, geo, persistent=True)
    _, src, _ = gen.generate()
    assert gen.tmem and gen.U == 6
    assert src.count("sf_tmem_alloc(") == 1 and src.count("sf_tmem_dealloc(") == 1
    assert src.index("sf_tmem_alloc(") < src.index("while (item <") < src.index("sf_tmem_dealloc(")
    # per unrolled step and field: one x8 + one x4 store and load of the 12 words; fast and boundary copies
    assert src.count("sf_tmem_st8(") == src.count("sf_tmem_ld8(") == 2 * 6 * 4
    assert src.count("sf_tmem_st4(") == src.count("sf_tmem_ld4(") == 2 * 6 * 4
    assert src.count("sf_tmem_wait_ld();") == 2 * 6 * 4
    # the switch off: the pass is what it was
    off = lower_stream.StreamKernelGen(prog, ops, ana, lower_stream.Geometry(ana, 4, 3, 24, 1, 5, 16),
                                       persistent=True).generate()[1]
    assert "sf_tmem" not in off


def _streamed(prog, **opts):
    from stencilflow_b200 import planner
    plan = planner.plan_program(prog, planner.PlanOptions(**opts) if opts else None)
    return [l for l in plan.lowered.launches if l.family == "streamed"]


def test_tmem_knob_reaches_the_generator():
    """diamond3d sits far below the register limit: tmem=1 keeps its planes in registers, tmem=2 parks them all the
    same, tmem=0 never parks; on the Jacobi-3D pass of config 1 (at its register limit) only tmem=0 keeps them."""
    geo = dict(max_depth=4, rows_per_thread=4, warps=8, threads_per_row=32, prefetch=2, sync="cta")
    prog = _program("diamond3d_12x10x16")
    assert [l.info["tmem"] for l in _streamed(prog, tmem=2, **geo)] == [{"a": 2, "r": 2}]
    assert [l.info["tmem_store"] for l in _streamed(prog, tmem=2, **geo)] == [{"a": 2, "r": -2}]
    assert [l.info["tmem"] for l in _streamed(prog, tmem=1, **geo)] == [{}]
    assert [l.info["tmem"] for l in _streamed(prog, tmem=0, **geo)] == [{}]
    # the register estimate, not the knob, decides at 1: 12 warps x 3 rows of config 1 parks, with the mbarriers
    config1 = dict(max_depth=4, rows_per_thread=3, warps=12, prefetch=5)
    prog = _program("ref_jacobi3d_32x32x32_8itr_8vec")
    on = _streamed(prog, tmem=1, **config1)
    assert [l.info["tmem"] for l in on] == [{"a": 2, "b0": 2, "b1": 2, "b2": 2}, {"b3": 2, "b4": 2, "b5": 2, "b6": 2}]
    assert all(l.info["sync"] == "flags" for l in on)
    assert not any(l.info["tmem"] for l in _streamed(prog, tmem=0, **config1))


def test_tmem_knob_from_the_environment(monkeypatch):
    from stencilflow_b200.planner import PlanOptions
    for value in ("0", "1", "2"):
        monkeypatch.setenv("SFB200_TMEM", value)
        assert PlanOptions().tmem == int(value) and not PlanOptions().is_default
    monkeypatch.delenv("SFB200_TMEM")
    assert PlanOptions().tmem == 1


@pytest.mark.parametrize("index,parked", [(1, True), (2, False), (3, False), (4, True)])
def test_default_plans_of_the_baseline_configs(monkeypatch, index, parked):
    """The cost model's policy: the Jacobi-3D passes of configs 1 and 4 park their planes and synchronise by
    per-field mbarriers; hdiff (config 2) and the 2-D chain (config 3) keep every plane in registers."""
    from stencilflow_b200 import programs
    from stencilflow_b200.planner import PlanOptions
    for knob in PlanOptions.KNOBS + ("SFB200_TUNED", "SFB200_PERSISTENT"):
        monkeypatch.delenv(knob, raising=False)
    name, prog, _ = programs.baseline_config(index)
    streamed = _streamed(_program_at(programs.write_program(prog, name)))
    assert streamed
    if parked:
        assert all(l.info["tmem"] and l.info["sync"] == "flags" for l in streamed)
    else:
        assert not any(l.info["tmem"] for l in streamed)


def test_gpu_matrix_covers_every_parking_shape(monkeypatch):
    """The GPU matrix of ``test_tmem_gpu.py``, lowered here: every entry parks what it says it parks, and together the
    entries reach every branch of the generator's parking code -- a slot parked at the start of the step (-2) and
    after an operator (>= 0), an age-3 slot, two fields parked at one point, float32 and float64, the chunk grid and
    persistent CTAs, and each synchronisation scheme.  Pruning the matrix must not drop one of them unnoticed."""
    import test_tmem_gpu as gm
    seen = set()
    for name, opts, env, slots in gm.MATRIX:
        for knob in ("SFB200_PERSISTENT", "SFB200_HALO_SKIP", "SFB200_SPLITLOOP"):
            monkeypatch.delenv(knob, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        prog = _program_at(gm.case_path(name))
        assert [l.info["tmem"] for l in _streamed(prog, tmem=0, **opts)] == [{}] * len(slots), (name, opts, env)
        on = _streamed(prog, tmem=2, **opts)
        assert [l.info["tmem"] for l in on] == slots, (name, opts, env)
        dtype = prog.ops[0].data_type.name
        for l in on:
            info = l.info
            if not info["tmem"]:
                continue
            points = list(info["tmem_store"].values())
            seen.update(("store", "start" if k == -2 else ("input" if k == -1 else "op")) for k in points)
            seen.update(("age", a) for a in info["tmem"].values())
            if len(points) > len(set(points)):
                seen.add("shared store point")
            seen.add(dtype)
            seen.add("persistent" if info["persistent"] else "chunk grid")
            seen.add(info["sync"])
            if info["direct"]:
                seen.add("direct")
            if info["halo_skip"][2] < len(l.ops):
                seen.add("halo warps")
    need = {("store", "start"), ("store", "op"), ("age", 1), ("age", 2), ("age", 3), "shared store point",
            "float32", "float64", "persistent", "chunk grid", "cta", "pair", "flags", "halves", "direct", "halo warps"}
    assert need <= seen, sorted(map(str, need - seen))


def test_chunk_grid_allocates_after_its_early_return(monkeypatch):
    """A CTA of the one-per-(tile, chunk) grid whose chunk is empty leaves before it allocates tensor memory; every
    other one frees its columns once, at the end."""
    from stencilflow_b200 import lower_stream
    monkeypatch.setenv("SFB200_PERSISTENT", "0")
    prog = _config1()
    ops = list(prog.ops)[:4]
    ana = _analysis(prog, ops)
    geo = lower_stream.Geometry(ana, 4, 3, 24, 1, 5, 16, "flags", tmem=True)
    gen = lower_stream.StreamKernelGen(prog, ops, ana, geo)
    _, src, _ = gen.generate()
    assert gen.tmem and not gen.persistent
    assert src.count("sf_tmem_alloc(") == 1 and src.count("sf_tmem_dealloc(") == 1
    assert src.index("if (c_begin >= c_end) return;") < src.index("sf_tmem_alloc(") < src.index("sf_tmem_dealloc(")
    assert "return;" not in src[src.index("sf_tmem_alloc("):]

"""Tensor-memory window slots of the fused 3-D pass (no GPU): which slots qualify, what the register estimate
and the shared-memory budget make of them, and what the generator emits."""
import pytest

from conftest import program_path


def _program(name):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    return make_program(KernelChainGraph(program_path(name)))


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

"""Host-side planning decisions (no GPU): the plans the BASELINE configs get, the options that reach
the generator, the chunking that fills every CTA slot of an SM."""
import os

import pytest

from conftest import program_path


def _program(index, variant=None):
    import bench
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    bench.VARIANT = variant
    try:
        name, prog, _ = bench.build_config(index)
    finally:
        bench.VARIANT = None
    return CudaProgram(programs.write_program(prog, name), allocate=False), prog


def test_config1_plan(native_lib):
    p, prog = _program(1)
    launches = p.lowered.launches
    assert [len(l.ops) for l in launches] == [4, 4] and all(l.family == "streamed" for l in launches)
    info = launches[0].info
    assert info["tile"] == [72, 64] and info["R"] == 3 and info["prefetch"] == 5 and info["unroll"] == 6
    assert launches[0].block == (384, 1, 1) and launches[0].smem <= 227 * 1024
    # persistent CTAs, one per SM, fetching items from a shared list: two waves of whole tiles, the 66
    # domain-edge tiles (slower: boundary code in every step) first, then the 8 tiles that do not fill a wave
    # in halving plane ranges so that the CTAs finish together
    assert info["persistent"] and info["tiles"] == 19 * 16
    assert launches[0].grid_fn(0, 1024) == (148, 1, 1)
    items = info["work_items_fn"](0, 1024)
    whole = items[:296]
    assert all((p0, p1) == (0, 1024) for _, p0, p1 in whole) and len({t for t, _, _ in whole}) == 296
    edge = {t for t in range(304) if t % 19 in (0, 18) or t // 19 in (0, 15)}
    assert {t for t, _, _ in whole[:len(edge)]} == edge
    rest = items[296:]
    assert len({t for t, _, _ in rest}) == 8 and not ({t for t, _, _ in rest} & {t for t, _, _ in whole})
    lengths = [p1 - p0 for _, p0, p1 in rest]
    assert lengths == sorted(lengths, reverse=True) and lengths[-1] <= 32
    for t in {t for t, _, _ in rest}:
        covered = sorted((p0, p1) for tt, p0, p1 in rest if tt == t)
        assert covered[0][0] == 0 and covered[-1][1] == 1024 and all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
    steps = sum(p1 - p0 + info["stream_overhead_planes"] for _, p0, p1 in items) / 148.0
    assert steps <= 1.02 * (19 * 16 * 1024 / 148.0)
    table = info["work_fn"](0, 1024)
    assert table[:3] == [0, 0, len(items)] and table[3:9] == [items[0][0], 0, 1024, items[1][0], 0, 1024]
    # algorithmic bytes of a pass: the field in, the field out
    assert launches[0].reads == ["a"] and launches[0].writes == ["b3"]


def test_config1_halving_list(native_lib, monkeypatch):
    """SFB200_SCHED=halving: the list the longest-first one replaced -- one wave of whole tiles (neighbours in
    lockstep), then the other 156 tiles in rounds of plane ranges that halve, 512, 256, ... 32."""
    monkeypatch.setenv("SFB200_SCHED", "halving")
    p, prog = _program(1)
    info = p.lowered.launches[0].info
    items = info["work_items_fn"](0, 1024)
    assert items[:148] == [(t, 0, 1024) for t in range(148)]
    rest = items[148:]
    assert {t for t, _, _ in rest} == set(range(148, 304))
    assert rest[:156] == [(t, 0, 512) for t in range(148, 304)]          # tile-minor: neighbours side by side
    lengths = [p1 - p0 for _, p0, p1 in rest]
    assert lengths == sorted(lengths, reverse=True) and lengths[-1] == 32
    for t in range(148, 304):
        covered = sorted((p0, p1) for tt, p0, p1 in rest if tt == t)
        assert covered[0][0] == 0 and covered[-1][1] == 1024 and all(a[1] == b[0] for a, b in zip(covered, covered[1:]))


@pytest.mark.parametrize("index", [1, 2, 3])
def test_cost_model_alone_finds_the_measured_plans(native_lib, monkeypatch, index):
    """SFB200_TUNED=0: without the table of measured plans the planner's cost model arrives at the same
    kernels for the three benchmark programs (the table is a record of measurements, not what the choice rests on)."""
    tuned = _program(index)[0]
    monkeypatch.setenv("SFB200_TUNED", "0")
    model = _program(index)[0]
    assert [l.kernel for l in model.lowered.launches] == [l.kernel for l in tuned.lowered.launches]
    assert [l.info["tile"] for l in model.lowered.launches] == [l.info["tile"] for l in tuned.lowered.launches]


def test_launch_bound_grids_are_not_fused(native_lib, tmp_path):
    """The latency terms of the cost model: on 32^3 ... 64^3 an 8-operator chain is eight one-operator launches
    (replayed through a CUDA graph), from 96^3 on it is fused passes (profiles/r02b_small_grid_sizes.txt)."""
    import json
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    for n, fused in ((32, False), (64, False), (96, True), (256, True)):
        path = tmp_path / "chain_{}.json".format(n)
        path.write_text(json.dumps(programs.jacobi3d_chain([n, n, n], 8)))
        p = CudaProgram(str(path), allocate=False)
        families = [l.family for l in p.lowered.launches]
        assert (families == ["streamed", "streamed"]) if fused else (families == ["general"] * 8), (n, families)


def test_pipelined_call_pieces_are_short_at_both_ends():
    """The overlapped host-array call: short pieces at both ends (what cannot overlap is the first upload and the
    last download), equal pieces in between, every plane exactly once."""
    from stencilflow_b200.cuda_program import CudaProgram
    for (n0, n1, pieces, reach) in [(0, 1024, 16, 4), (0, 32768, 16, 8), (100, 612, 8, 2), (0, 80, 16, 1), (0, 2048, 32, 4)]:
        ends = CudaProgram._piece_ends(n0, n1, pieces, reach)
        sizes = [b - a for a, b in zip([n0] + ends[:-1], ends)]
        assert ends[-1] == n1 and all(s_ > 0 for s_ in sizes) and ends == sorted(ends)
        if (n1 - n0) // pieces > 8 * reach:
            assert sizes[0] == max(4 * reach, 8) == sizes[-1] and sizes[0] < max(sizes)
            assert sizes[1] == 2 * sizes[0] == sizes[-2] and sizes == sizes[::-1][:len(sizes)] or sum(sizes) == n1 - n0
            assert sum(1 for s_ in sizes if s_ >= max(sizes) - 1) >= pieces // 2
    os.environ["SFB200_PIPELINE_RAMP"] = "0"
    try:
        assert CudaProgram._piece_ends(0, 1024, 16, 4) == [64 * (s_ + 1) for s_ in range(16)]
    finally:
        del os.environ["SFB200_PIPELINE_RAMP"]


def test_config3_plan_uses_small_independent_ctas(native_lib, monkeypatch):
    p, prog = _program(3)
    launches = p.lowered.launches
    assert [len(l.ops) for l in launches] == [8, 8]
    l = launches[0]
    # one-warp CTAs, eight of them per SM (255 registers each), each with its own TMA ring and barrier
    assert l.block == (32, 1, 1) and l.info["tile"] == [1, 128] and l.info["prefetch"] == 5
    # 293 column tiles on 8 x 148 CTA slots: fewer tiles than slots, so the plain (tile, chunk) grid is used
    assert not l.info["persistent"] and l.info["tiles"] == 293
    gx, gy, gz = l.grid_fn(0, 32768)
    assert gx == 293 and gy == 1
    # many short chunks (at most 32 x the 16 warm-up rows each: measured 4.7 % faster than the few long chunks
    # that minimise waves x (rows + warm-up)), the last wave of CTAs nearly full
    waves = gx * gz / (8 * 148.0)
    assert waves >= 12 and (waves - int(waves) > 0.8 or waves == int(waves))
    assert l.info["chunk_fn"](0, 32768) <= 32 * l.info["stream_overhead_planes"]
    assert l.info["stream_overhead_planes"] * gz <= 0.04 * 32768
    # ... unless persistent CTAs are forced: every tile cut into row ranges, long ones first
    monkeypatch.setenv("SFB200_PERSISTENT", "1")
    p, prog = _program(3)
    l = p.lowered.launches[0]
    items = l.info["work_items_fn"](0, 32768, 8 * 148)
    assert l.info["persistent"] and l.grid_fn(0, 32768, 8 * 148) == (min(8 * 148, len(items)), 1, 1)
    assert [t for t, _, _ in items[:293]] == list(range(293))          # tile-minor: neighbours side by side
    rows = sorted((p0, p1) for (t, p0, p1) in items if t == 5)
    assert rows[0][0] == 0 and rows[-1][1] == 32768 and all(a[1] == b[0] for a, b in zip(rows, rows[1:]))
    overhead = l.info["stream_overhead_planes"]
    assert min(p1 - p0 for p0, p1 in rows) >= 4 * overhead


def test_one_cta_per_tile_chunk_grid_still_available(native_lib, monkeypatch):
    monkeypatch.setenv("SFB200_PERSISTENT", "0")
    p, prog = _program(1)
    l = p.lowered.launches[0]
    assert not l.info["persistent"] and ("chunk",) in l.args
    gx, gy, gz = l.grid_fn(0, 1024)
    assert (gx, gy) == (19, 16) and gx * gy * gz >= 4 * 148


@pytest.mark.parametrize("sched", ["lpt", "rows", "halving"])
def test_schedule_work_covers_every_plane_once(monkeypatch, sched):
    from stencilflow_b200.lower_stream import schedule_work, pack_work_table
    monkeypatch.setenv("SFB200_SCHED", sched)
    for (tiles, planes, slots, ov) in [(304, 1024, 148, 8), (1184, 256, 148, 8), (150, 1024, 148, 8), (1, 32, 148, 8),
                                       (24, 1024, 148, 5), (137, 32768, 592, 16), (3, 7, 148, 2), (600, 64, 148, 8),
                                       (304, 64, 148, 8), (2, 1024, 148, 8), (1184, 2048, 148, 8), (296, 1024, 148, 8),
                                       (297, 40, 148, 8)]:
        # (domain-edge tiles as the lowering passes them: a frame around a 19-wide grid of tiles)
        edge = {t for t in range(tiles) if t % 19 in (0, 18) or t < 19 or t >= tiles - 19}
        items = schedule_work(tiles, planes, slots, ov, edge_tiles=edge)
        seen = {}
        for (t, p0, p1) in items:
            assert 0 <= t < tiles and 0 <= p0 < p1 <= planes
            seen.setdefault(t, []).append((p0, p1))
        assert sorted(seen) == list(range(tiles))
        for t, ranges in seen.items():
            ranges.sort()
            assert ranges[0][0] == 0 and ranges[-1][1] == planes
            assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        # longest items first: what is fetched late is short
        lengths = [p1 - p0 for _, p0, p1 in items]
        assert lengths[0] == max(lengths)
        # the warm-up planes every item re-streams stay a small part of a big pass
        if tiles * planes >= 64 * slots * ov:
            assert sum(p1 - p0 + ov for _, p0, p1 in items) <= 1.06 * tiles * planes
        table = pack_work_table(items)
        assert table[:3] == [0, 0, len(items)] and len(table) == 3 + 3 * len(items)
    # exactly 8 tiles per SM (config 4 on 8 GPUs): whole tiles only, nothing is cut
    assert schedule_work(1184, 256, 148, 8) == [(t, 0, 256) for t in range(1184)]
    # a tiny grid is cut as finely as its single tile allows: launch latency, not warm-up, is what counts
    assert len(schedule_work(1, 32, 148, 8)) == 32


def test_cost_model_picks_small_ctas_and_depth_for_untuned_2d(native_lib):
    p, prog = _program(3, "w1d")                      # not in the table of measured plans
    launches = p.lowered.launches
    assert [len(l.ops) for l in launches] == [8, 8]
    assert launches[0].block == (32, 1, 1) and launches[0].info["prefetch"] == 5     # one-warp CTAs, eight per SM
    assert "w" in launches[0].reads                   # the 1-D weight is read by the fused pass itself


def test_direct_rows_option_reaches_the_generator(native_lib):
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    path = program_path("ref_jacobi3d_32x32x32_8itr_8vec")
    on = CudaProgram(path, allocate=False, plan_options=PlanOptions(max_depth=4, rows_per_thread=4, warps=8,
                                                                     threads_per_row=32, prefetch=4, direct=1))
    off = CudaProgram(path, allocate=False, plan_options=PlanOptions(max_depth=4, rows_per_thread=4, warps=8,
                                                                      threads_per_row=32, prefetch=4))
    assert on.lowered.launches[0].info["direct"] == ["a"] and off.lowered.launches[0].info["direct"] == []
    # no exchange ring for the input, one more TMA slot instead
    src_on = on.lowered.kernels[on.lowered.launches[0].kernel].source
    src_off = off.lowered.kernels[off.lowered.launches[0].kernel].source
    assert "xrow_f0" not in src_on and "xrow_f0" in src_off
    # a non-zero boundary value needs the fix-up in registers: the option leaves that input on the ring
    keep = CudaProgram(program_path("jacobi3d_16x24x32_5itr_const1"), allocate=False,
                       plan_options=PlanOptions(max_depth=4, rows_per_thread=4, warps=8, threads_per_row=32,
                                                prefetch=4, direct=1))
    assert keep.lowered.launches[0].info["direct"] == []


def test_environment_knobs(monkeypatch):
    from stencilflow_b200.planner import PlanOptions
    for k in PlanOptions.KNOBS:
        monkeypatch.delenv(k, raising=False)
    assert PlanOptions().is_default
    monkeypatch.setenv("SFB200_DIRECT", "1")
    monkeypatch.setenv("SFB200_SYNC", "pair")
    o = PlanOptions()
    assert o.direct == 1 and o.sync == "pair" and not o.is_default
    assert PlanOptions(direct=0).direct == 0


def test_reference_arm_line(monkeypatch):
    """`bench.py --impl reference`: one JSON line with the contract's keys, timed on all host threads
    even when the launcher exports OMP_NUM_THREADS=1 (torchrun does), the thread count taken from the
    OpenMP runtime itself."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    env = dict(os.environ, OMP_NUM_THREADS="1")
    env.pop("SFB200_REF_THREADS", None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "0",
                          "--steps", "3", "--warmup", "1"], stdout=subprocess.PIPE, text=True, env=env, timeout=300,
                         check=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "stencil_cell_updates_per_s"
    assert line["unit"] == "cell-updates/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["ms_per_step"] > 0 and "32x32x32" in line["config"]["workload"]
    # exactly the requested number of timed executions; the same config keys as the GPU arm prints
    assert line["steps"] == 3 and line["warmup"] == 1
    assert set(line["config"]) == {"workload", "per_gpu", "l2", "input"}


def test_bench_dump_outputs_writes_a_fixed_sample(tmp_path):
    """``bench.py --dump-outputs``: a small output is written whole, a large one as the same seeded sample
    on every run, all files within the size budget; the undefined -halo border is left out."""
    import types
    import numpy as np
    import bench
    fields = {"small": np.arange(6 * 7 * 8, dtype=np.float64).reshape(6, 7, 8),
              "large": np.full((68, 512, 260), np.nan, np.float32)}
    fields["large"][2:-2, 2:-2, 2:-2] = np.random.default_rng(0).random((64, 508, 256), np.float32)
    fake = types.SimpleNamespace(program=types.SimpleNamespace(outputs=list(fields)),
                                 download=lambda name: fields[name].copy())
    for run in ("a", "b"):
        bench.dump_outputs(fake, str(tmp_path / run), halo=2)
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), fields["small"][2:-2, 2:-2, 2:-2])
    large = np.load(tmp_path / "a" / "large.npy")
    assert large.dtype == np.float32 and large.ndim == 1 and large.size > 1000000
    assert not np.isnan(large).any()
    assert np.array_equal(large, np.load(tmp_path / "b" / "large.npy"))
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 << 20


def test_choose_chunk_balances_waves_and_warmup():
    from stencilflow_b200.lower_stream import choose_chunk
    # 304 tiles of config 1, 8 warm-up planes per chunk, one CTA per SM
    ci = choose_chunk(1024, 304, 8, sms=148)

    def cost(c):                                  # rounds of CTAs x planes each CTA streams
        return -(-(304 * -(-1024 // c)) // 148) * (c + 8)
    assert cost(ci) == min(cost(-(-1024 // n)) for n in range(1, 65)) and 8.0 / ci < 0.08
    # a single tile column must be cut into many chunks to occupy the machine at all
    ci = choose_chunk(32768, 1, 16, sms=148)
    assert -(-32768 // ci) >= 60
    # more resident CTAs per SM -> more, shorter chunks
    assert choose_chunk(32768, 137, 16, sms=4 * 148) < choose_chunk(32768, 137, 16, sms=148)


@pytest.mark.parametrize("name,depth,expect", [
    ("ref_jacobi3d_32x32x32_8itr_8vec", 4, (4, 8)),      # two passes of four: 4 per pass, 8 in total
    ("ref_jacobi3d_32x32x32_8itr_8vec", 2, (2, 8)),
    ("ref_jacobi3d_32x32x32_8itr_8vec", 8, (8, 8)),
    ("hdiff_24x28x16", 4, (2, 2)),                        # lap -> flx/fly -> out reaches 2 planes along i
])
def test_halo_depth_and_total_reach(native_lib, name, depth, expect):
    from stencilflow_b200 import distributed
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    p = CudaProgram(program_path(name), allocate=False, plan_options=PlanOptions(max_depth=depth))
    assert (distributed.halo_depth(p.lowered), distributed.total_reach(p.lowered)) == expect


def test_halo_schedule_of_a_two_pass_chain(native_lib):
    from stencilflow_b200 import distributed
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    p = CudaProgram(program_path("ref_jacobi3d_32x32x32_8itr_8vec"), allocate=False,
                    plan_options=PlanOptions(max_depth=4))
    middle = distributed.Slab(1, 4, 32, 4)
    sends = distributed.halo_schedule(p.lowered, middle)
    # only the first pass's result crosses slab boundaries: 4 planes up, 4 planes down
    assert sorted((s.launch, s.field, s.peer, s.src_end - s.src_begin) for s in sends) == \
        [(0, "b3", 0, 4), (0, "b3", 2, 4)]
    assert distributed.halo_schedule(p.lowered, distributed.Slab(0, 1, 32, 4)) == []


def test_partition_cache_distinguishes_source_type(native_lib, tmp_path):
    """Two chains with identical taps but sources of different type: float32 operators on a float32
    field stream, the same operators on a float64 field cannot (mixed types) -- the cost cache of the
    partition must not carry the first answer over to the second (either order)."""
    import json
    from stencilflow_b200.cuda_program import CudaProgram

    def chain(src, names):
        out, prev = {}, src
        for n in names:
            out[n] = {"data_type": "float32", "boundary_conditions": {prev: {"type": "constant", "value": 0.0}},
                      "computation_string": "{n} = 0.25 * ({p}[i,j,k-1] + {p}[i,j,k+1] + {p}[i-1,j,k] + {p}[i,j+1,k])".format(n=n, p=prev)}
            prev = n
        return out

    for order in ((("a", "float32"), ("b", "float64")), (("b", "float64"), ("a", "float32"))):
        prog = {"dimensions": [96, 128, 256], "outputs": [], "inputs": {}, "program": {}}
        for k, (src, dt) in enumerate(order):
            prog["inputs"][src] = {"data": "constant:1.0", "data_type": dt}
            names = ["o{}_{}".format(src, s) for s in range(3)]
            prog["program"].update(chain(src, names))
            prog["outputs"].append(names[-1])
        path = tmp_path / "mixed_{}.json".format(order[0][0])
        path.write_text(json.dumps(prog))
        p = CudaProgram(str(path), allocate=False)            # must plan without raising in either order
        fam = {op: l.family for l in p.lowered.launches for op in l.ops}
        group = {op: tuple(l.ops) for l in p.lowered.launches for op in l.ops}
        # the float32 chain on the float32 field streams (its first stage may be cheaper as a one-operator
        # launch on a grid this small: a streamed kernel costs a few microseconds before its first plane) ...
        assert all(fam["oa_{}".format(k)] == "streamed" for k in (1, 2)), (fam, group)
        # ... the operator reading the float64 field into a float32 result cannot (mixed types)
        assert fam["ob_0"] == "general", (fam, group)

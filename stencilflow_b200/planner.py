"""Fusion-depth and tile planner: decides how the operator DAG is cut into passes over HBM.

This replaces the reference's buffer-placement optimizer (``stencilflow/optimizer.py:73-307``), which
greedily moves FPGA delay/window buffers between fast (on-chip) and slow (off-chip) memory under a
size or communication-volume bound.  On a GPU the same trade-off reads: a field that stays *inside* a
pass lives in registers/shared memory (fast memory) and costs no HBM traffic; a field that crosses a
pass boundary is written to and re-read from HBM (slow memory).  The planner therefore

1. walks the operators in topological order and grows a *pass* (fusion group) while the group is
   streamable (see :mod:`lower_stream` for the conditions), its fusion depth stays within
   ``max_depth`` and its tile fits the shared-memory/register budget (227 KB per CTA, 64 K registers
   per SM);
2. lowers each pass with the streamed template, or -- for operators the template cannot express
   (copy boundaries, far taps, lower-dimensional array inputs, mixed boundary values ...) -- with the
   general one-operator kernel;
3. assigns HBM storage to the fields that cross pass boundaries, reusing the storage of dead
   intermediates (the reference keeps every transient alive, ``stencilflow/sdfg_generator.py:626-630``;
   results are identical, the footprint is what makes 2048^3 x 64 operators fit).

``Plan.describe()`` is the inspectable record of these decisions (written to ``plan.json`` next to
the generated source).
"""

import hashlib
import json
import os
from typing import Dict, List, Optional

from . import lower_cuda
from .stencil_op import StencilProgram


# default of PlanOptions.tmem (SFB200_TMEM): park window planes in tensor memory where a 3-D pass needs the registers
TMEM_DEFAULT = "1"
TUNED_PLANS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tuned_plans.json")


def structure_key(program: StencilProgram) -> str:
    """Hash of the operator structure that determines the best plan, independent of names, extents
    and chain length: the *set* of distinct operator signatures, an operator's signature being its
    type, its boundary handling and its taps with each source named relative to the operator (the
    n-th operator before it, or the n-th program input).  An 8- and a 64-stage chain of the same
    stencil share a key; ``lookup_tuned`` then picks the entry with the closest extents."""
    op_index = {op.name: n for n, op in enumerate(program.ops)}
    inputs = [name for name, f in program.fields.items() if f.kind == "input"]

    def rel(field, k):
        if field in op_index:
            return "op-{}".format(k - op_index[field])
        return "in{}".format(inputs.index(field)) if field in inputs else field

    sigs = set()
    for k, op in enumerate(program.ops):
        taps = sorted((rel(f, k), tuple(map(tuple, op.offsets3(f)))) for f in op.accesses)
        bcs = sorted((rel(f, k), bc.get("btype"), repr(bc.get("value")))
                     for f, bc in op.boundary_conditions.items() if f in op.accesses)
        sigs.add(json.dumps([op.data_type.name, taps, bcs, len(op.statements)], default=str))
    text = json.dumps([len(program.shape), sorted(sigs)])
    return hashlib.sha1(text.encode()).hexdigest()[:16]


def lookup_tuned(program: StencilProgram, table=None):
    """Entry of the measured-plan table for ``program``: same operator structure, and the extents
    closest (in log distance) among the entries whose innermost dimension is in the same class
    (narrow / wide) and whose cell count is within 64x.  None if there is none."""
    import math
    table = load_tuned() if table is None else table
    entries = table.get(structure_key(program))
    if not entries:
        return None
    shape = list(program.shape)
    best = None
    for entry in entries:
        other = entry.get("shape")
        if not other or len(other) != len(shape) or (other[-1] < 128) != (shape[-1] < 128):
            continue
        dist = sum(abs(math.log2(a / float(b))) for a, b in zip(shape, other))
        if dist > 6.0:
            continue
        if best is None or dist < best[0]:
            best = (dist, entry)
    return best[1] if best else None


def load_tuned():
    """The table ``scripts/tune.py`` measures on a B200: structure key -> plan options."""
    try:
        with open(TUNED_PLANS) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


class PlanOptions:
    """Knobs, all overridable through ``SFB200_*`` environment variables.  When neither the caller
    nor the environment sets any of them, ``plan_program`` looks the program up in the table of
    measured plans (``tuned_plans.json``) before falling back on the cost model."""

    KNOBS = ("SFB200_FUSE", "SFB200_MAX_DEPTH", "SFB200_ROWS", "SFB200_WARPS", "SFB200_CHUNK", "SFB200_PREFETCH",
             "SFB200_VEC", "SFB200_KS", "SFB200_SYNC", "SFB200_DIRECT",
             "SFB200_TMEM")

    def __init__(self, fuse=None, max_depth=None, rows_per_thread=None, warps=None, chunk=None,
                 prefetch=None, vector=None, threads_per_row=None, sync=None, direct=None, tmem=None,
                 peer_push=None, cluster=None, unaligned=None):
        env = os.environ
        self.is_default = (all(v is None for v in (fuse, max_depth, rows_per_thread, warps, chunk, prefetch, vector,
                                                   threads_per_row, sync, direct, tmem))
                           and not any(k in env for k in self.KNOBS) and env.get("SFB200_TUNED", "1") != "0")
        self.vector = int(env.get("SFB200_VEC", "0")) if vector is None else vector
        self.threads_per_row = int(env.get("SFB200_KS", "0")) if threads_per_row is None else threads_per_row
        self.fuse = (env.get("SFB200_FUSE", "1") != "0") if fuse is None else fuse
        self.max_depth = int(env.get("SFB200_MAX_DEPTH", "0")) if max_depth is None else max_depth
        self.rows_per_thread = int(env.get("SFB200_ROWS", "0")) if rows_per_thread is None else rows_per_thread
        self.warps = int(env.get("SFB200_WARPS", "0")) if warps is None else warps
        self.chunk = int(env.get("SFB200_CHUNK", "0")) if chunk is None else chunk
        self.prefetch = int(env.get("SFB200_PREFETCH", "0")) if prefetch is None else prefetch
        self.sync = env.get("SFB200_SYNC", "") if sync is None else sync
        # 1: neighbour rows of a streamed *input* field are read straight from its TMA ring (which then
        # keeps a plane one step longer) instead of being re-published through an exchange ring
        self.direct = int(env.get("SFB200_DIRECT", "0")) if direct is None else int(direct)
        # 1: 3-D passes with one CTA per SM that sit at their register limit park the oldest plane of a window in
        # tensor memory between its last use as a centre plane and its use as an own-cell operand; 2: park every
        # slot that qualifies, whatever the register estimate (tests); 0: never
        self.tmem = int(env.get("SFB200_TMEM", TMEM_DEFAULT)) if tmem is None else int(tmem)
        # 1: a program whose fields fit the distributed shared memory of one 8-CTA cluster runs as one launch of
        # the cluster family (lower_cluster); 0: never.  Like ``peer_push`` not a tuning knob: it does not take
        # part in ``is_default`` and survives the replacement of the options by a measured plan.  Ignored with
        # fuse=False and in slab mode.
        self.cluster = int(env.get("SFB200_CLUSTER", "0")) if cluster is None else int(cluster)
        # 1: groups whose innermost row is not a multiple of 16 bytes stream too: the threads copy their input cells
        # into the shared-memory ring with cp.async (a tiled TMA map needs 16-byte row strides), and results leave by
        # single-cell stores (lower_stream).  0: such groups run as one-operator kernels.  Programs with aligned rows
        # get the same kernels either way.  Like ``cluster`` not a tuning knob; ignored with fuse=False and in slab mode.
        self.unaligned = int(env.get("SFB200_UNALIGNED", "0")) if unaligned is None else int(unaligned)
        # slab mode (set by distributed.SlabProgram): streamed kernels store the edge planes of their
        # results straight into the neighbouring GPUs' halo planes.  Not a tuning knob: it does not
        # take part in ``is_default`` and survives the replacement of the options by a measured plan.
        self.peer_push = bool(peer_push)

    def as_dict(self):
        return {k: v for k, v in self.__dict__.items() if k != "is_default"}


def share_storage(steps, nbytes, own=()) -> Dict[str, int]:
    """field -> storage id for the fields written by ``steps``, a sequence of (reads, writes) in execution
    order.  The fields in ``own`` come first, each with storage of its own.  Every other field takes the
    storage of a field of the same byte size that no step at or after its own writer reads, else new
    storage."""
    last_read = {}
    for idx, (reads, writes) in enumerate(steps):
        for f in reads:
            last_read[f] = idx
    assign, next_id = {}, 0
    free_pool = []            # (nbytes, storage id)
    busy = []                 # (last read index, nbytes, storage id)
    for name in own:
        assign[name] = next_id
        next_id += 1
    for idx, (reads, writes) in enumerate(steps):
        still = []
        for (lr, nb, sid) in busy:
            if lr < idx:
                free_pool.append((nb, sid))
            else:
                still.append((lr, nb, sid))
        busy = still
        for f in writes:
            if f in assign:
                continue
            nb = nbytes[f]
            sid = None
            for k, (pnb, psid) in enumerate(free_pool):
                if pnb == nb:
                    sid = psid
                    free_pool.pop(k)
                    break
            if sid is None:
                sid = next_id
                next_id += 1
            assign[f] = sid
            busy.append((last_read.get(f, idx), nb, sid))
    return assign


class Plan:
    def __init__(self, program: StencilProgram, lowered, passes, options):
        self.program = program
        self.lowered = lowered
        self.passes = passes          # list of dicts: {"ops": [...], "family": ..., ...}
        self.options = options

    def materialized_fields(self) -> List[str]:
        names = []
        for l in self.lowered.launches:
            for f in list(l.reads) + list(l.writes):
                if f not in names and not self.program.fields[f].is_scalar:
                    names.append(f)
        for name, f in self.program.fields.items():
            if f.kind in ("input", "output") and not f.is_scalar and name not in names:
                names.append(name)
        return names

    def buffer_assignment(self) -> Dict[str, int]:
        """field -> storage id.  Inputs and outputs own their storage; intermediates that cross
        pass boundaries share storage once dead (equal byte size only)."""
        fields = self.program.fields
        own = [name for name in self.materialized_fields() if fields[name].kind != "intermediate"]
        return share_storage([(l.reads, l.writes) for l in self.lowered.launches],
                             {name: f.nbytes for name, f in fields.items()}, own)

    def algorithmic_bytes(self) -> int:
        return self.lowered.algorithmic_bytes()

    def cell_updates(self) -> int:
        return len(self.program.ops) * self.program.cells

    def describe(self):
        fields = self.program.fields
        return {
            "program": self.program.name,
            "shape": list(self.program.shape),
            "operators": len(self.program.ops),
            "cell_updates": self.cell_updates(),
            "options": self.options.as_dict(),
            "tuned_from": getattr(self, "tuned_from", None),
            "passes": [
                {
                    "family": l.family, "kernel": l.kernel, "ops": l.ops, "reads": l.reads,
                    "writes": l.writes, "block": list(l.block), "smem": l.smem,
                    "algorithmic_bytes": sum(fields[f].nbytes for f in l.reads) +
                    sum(fields[f].nbytes for f in l.writes),
                    "info": {k: v for k, v in l.info.items() if not callable(v)},
                } for l in self.lowered.launches
            ],
            "algorithmic_bytes": self.algorithmic_bytes(),
            "storage": self.buffer_assignment(),
        }


def plan_program(program: StencilProgram, options: Optional[PlanOptions] = None,
                 specialize=None) -> Plan:
    options = options or PlanOptions()
    tuned_from = None
    if options.is_default:
        entry = lookup_tuned(program)
        if entry:
            options = PlanOptions(**dict(entry["options"], peer_push=options.peer_push, cluster=options.cluster,
                                         unaligned=options.unaligned))
            tuned_from = entry.get("measured")
    lowered = lower_cuda.LoweredProgram(program)
    passes = []
    groups = None
    if options.cluster and options.fuse and not options.peer_push:
        from . import lower_cluster
        layout = lower_cluster.ClusterLayout(program)
        if layout.fits:
            lower_cluster.lower_program_cluster(lowered, layout, specialize)
            plan = Plan(program, lowered, [{"family": "cluster", "ops": [op.name for op in program.ops]}], options)
            plan.tuned_from = tuned_from
            return plan
    if options.fuse:
        try:
            from . import lower_stream
        except ImportError:
            lower_stream = None
        if lower_stream is not None:
            groups = lower_stream.partition(program, options)
    if groups is None:
        groups = [("general", [op]) for op in program.ops]
    for family, ops in groups:
        if family == "general":
            for op in ops:
                lower_cuda.lower_general_op(lowered, op, specialize)
                passes.append({"family": "general", "ops": [op.name]})
        else:
            from . import lower_stream
            try:
                lower_stream.lower_group(lowered, ops, options, specialize)
                passes.append({"family": "streamed", "ops": [op.name for op in ops]})
            except lower_stream.NotStreamable:
                # the partition's estimate was wrong about this group: one-operator kernels always work
                for op in ops:
                    lower_cuda.lower_general_op(lowered, op, specialize)
                    passes.append({"family": "general", "ops": [op.name]})
    plan = Plan(program, lowered, passes, options)
    plan.tuned_from = tuned_from
    return plan

"""The ``cluster`` kernel family: a whole small program in one launch of one thread-block cluster.

Grids of a few thousand cells are bound by launch latency, not by any pipe (DESIGN §3.4).  When every
field the program keeps fits the distributed shared memory of one cluster of C <= 8 CTAs (the portable
cluster size), all operators run in one kernel:

* **Ownership.** The outermost dimension (i in 3-D, j in 2-D, k in 1-D) is cut into C contiguous
  ranges of P planes (rows, or k-cells that are a multiple of the widest vector), one per CTA.  A CTA
  holds its range of every field that lives in shared memory, at the same offset in every CTA.
* **Shared memory.** Full-dimensional inputs are copied from HBM into the owner's shared memory once, at
  kernel start.  Results read by a later operator stay in shared memory; slots are reused once a field is
  dead (:func:`planner.share_storage`).  Lower-dimensional and 0-D inputs are read as ``sf_general``
  reads them: global memory and kernel arguments.
* **Operators** run in topological order, each CTA computing its own cells, V consecutive k-cells per
  thread.  The per-cell code is :meth:`GeneralKernelGen.emit_cell` -- the same tap grouping, boundary
  selects, compute type, literals and statements -- so the results are bit-identical to the one-operator
  kernels.  Only the row source differs: a row of another CTA is addressed through ``mapa`` (distributed
  shared memory), a row of the thread's own range is a local shared-memory address.
* **Synchronisation.** A cluster barrier (release/acquire) goes before an operator that reads a field
  written, or writes a slot read or written, since the previous barrier; one more precedes the exit so
  that no CTA leaves while a peer still reads its shared memory.

The cluster size is compile-time (``__cluster_dims__``), so the launch is a plain ``cuLaunchKernel`` of
grid (C, 1, 1).
"""

import hashlib

from .lower_cuda import GeneralKernelGen, KernelSpec, LaunchSpec, ctype_of, vector_width

CLUSTER_MAX = 8                  # portable cluster size
SMEM_LIMIT = 227 * 1024          # dynamic shared memory a CTA may opt into on sm_100a
MAX_THREADS = 1024
MAX_ITEMS_PER_THREAD = 8         # V-cell items a thread computes per operator (48^3 Jacobi-3D: 3.4)
SLOT_ALIGN = 16

CLUSTER_PRELUDE = r"""
// ---- thread-block cluster / distributed shared memory (sm_90+) ----
__device__ __forceinline__ u32 sf_cluster_rank() {
    u32 r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// generic address of the same shared-memory variable in CTA `rank` of the cluster
template <typename T>
__device__ __forceinline__ const T* sf_cl_map(const T* p, u32 rank) {
    u64 r;
    asm("mapa.u64 %0, %1, %2;" : "=l"(r) : "l"(p), "r"(rank));
    return reinterpret_cast<const T*>(r);
}
// element k of a 1-D field cut into chunks of P cells, one per CTA (an out-of-range k is never dereferenced;
// it is clamped so that the address handed to mapa stays inside a slot)
template <typename T, int P, int C>
__device__ __forceinline__ const T* sf_cl_at(const T* slot, int k) {
    const int kc = min(max(k, 0), C * P - 1);
    const int o = kc / P;
    return sf_cl_map(slot + (kc - o * P), (u32)o);
}
// a 0-D input as the loop body sees it: opaque, so that nothing computed from it alone is hoisted out of the
// loop over a thread's cells (a product of two scalars computed once before the loop is rounded on its own,
// where the one-operator kernel contracts it into an FMA with the sum it belongs to)
__device__ __forceinline__ float sf_keep(float x) { asm volatile("" : "+f"(x)); return x; }
__device__ __forceinline__ double sf_keep(double x) { asm volatile("" : "+d"(x)); return x; }
__device__ __forceinline__ int sf_keep(int x) { asm volatile("" : "+r"(x)); return x; }
__device__ __forceinline__ unsigned sf_keep(unsigned x) { asm volatile("" : "+r"(x)); return x; }
__device__ __forceinline__ long long sf_keep(long long x) { asm volatile("" : "+l"(x)); return x; }
__device__ __forceinline__ unsigned long long sf_keep(unsigned long long x) { asm volatile("" : "+l"(x)); return x; }
template <typename T>
__device__ __forceinline__ T sf_keep(T x) { return (T)sf_keep((int)x); }
__device__ __forceinline__ void sf_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
"""


def _ceil(a, b):
    return -(-a // b)


class ClusterLayout:
    """Host-side plan of a cluster kernel: ownership, shared-memory slots, barriers and block size.
    ``fits`` is the capacity rule (checked before any code is generated)."""

    def __init__(self, program):
        from .planner import share_storage
        self.program = program
        fields = program.fields
        ops = program.ops
        self.outer = program.iterators[0]
        self.n = program.shape[0]
        self.vecs = [vector_width(program, op) for op in ops]
        unit = max(self.vecs) if len(program.shape) == 1 else 1
        units = self.n // unit
        c = min(CLUSTER_MAX, units)
        p_units = _ceil(units, c)
        self.C = _ceil(units, p_units)                   # fewer CTAs if the last ranges would be empty
        self.P = p_units * unit                          # planes / rows / k-cells per CTA
        self.plane = program.cells // self.n             # elements per index of the outermost dimension
        self.ranges = [[c * self.P, min(self.n, (c + 1) * self.P)] for c in range(self.C)]
        full = list(program.iterators)
        read_later = {f for op in ops for f in op.accesses}
        self.inputs = [name for name, f in fields.items()
                       if f.kind == "input" and not f.is_scalar and name in read_later]
        self.loaded = [name for name in self.inputs if fields[name].dims == full]
        self.smem = self.loaded + [op.name for op in ops if op.name in read_later]
        slot_bytes = {f: _ceil(self.P * self.plane * fields[f].data_type.bytes, SLOT_ALIGN) * SLOT_ALIGN
                      for f in self.smem}
        steps = [([], list(self.loaded))]
        steps += [([f for f in op.accesses if f in slot_bytes], [op.name] if op.name in slot_bytes else [])
                  for op in ops]
        sid = share_storage(steps, slot_bytes)
        offsets, total = {}, 0
        for s in sorted(set(sid.values())):
            offsets[s] = total
            total += next(slot_bytes[f] for f in sid if sid[f] == s)
        self.slot = {f: sid[f] for f in self.smem}
        self.offset = {f: offsets[sid[f]] for f in self.smem}
        self.smem_bytes = total
        # barriers: before op m when it reads a field written, or writes a slot read or written, since the last one
        self.barriers = []
        written, touched = set(self.loaded), set()
        for m, op in enumerate(ops):
            reads = [f for f in op.accesses if f in self.slot]
            mine = self.slot.get(op.name)
            if any(f in written for f in reads) or (mine is not None and (
                    mine in touched or mine in {self.slot[f] for f in written})):
                self.barriers.append(m)
                written, touched = set(), set()
            touched |= {self.slot[f] for f in reads}
            if mine is not None:
                written.add(op.name)
        items = max(_ceil(self.P * self.plane, v) for v in self.vecs)
        self.threads = min(MAX_THREADS, _ceil(items, 32) * 32)
        # capacity: the CTA's slots fit its shared memory, and its cells fit a few items per thread (a program that
        # keeps nothing in shared memory must not run a large grid on C SMs)
        self.fits = self.smem_bytes <= SMEM_LIMIT and items <= MAX_ITEMS_PER_THREAD * MAX_THREADS

    def describe(self):
        return {"cluster": self.C, "outer": self.outer, "planes_per_cta": self.P, "ranges": self.ranges,
                "slots": {f: [self.offset[f], self.slot[f]] for f in self.smem}, "barriers_before": self.barriers,
                "threads": self.threads}


class ClusterOpGen(GeneralKernelGen):
    """One operator's per-cell code inside the cluster kernel: rows of fields in shared memory come
    from the owning CTA; everything else is the general kernel's."""

    def __init__(self, op, program, layout, specialize=None):
        super().__init__(op, program, specialize)
        self.layout = layout
        self.slab_axis = None           # one cluster computes the whole domain

    def _row_pointer(self, field, di, dj, rid, base):
        lay = self.layout
        if field not in lay.slot:
            return super()._row_pointer(field, di, dj, rid, base)
        ft = ctype_of(self.program.fields[field].data_type)
        slot = "sm{}".format(lay.smem.index(field))
        NI, NJ, NK = self.n3
        if lay.outer == "k":
            return "  const {}* __restrict__ p{} = {};".format(ft, rid, slot)
        if lay.outer == "i":
            pos, off, rest = "i", di, " + (j + ({})) * {}".format(dj, NK)
        else:
            pos, off, rest = "j", dj, ""
        if not off:
            return "  const {}* __restrict__ p{} = {} + ({} - lo) * {}{};".format(ft, rid, slot, pos, lay.plane, rest)
        # a masked row is never read, but the address handed to mapa stays inside the owner's slot: the row
        # falls back to the thread's own (i, j)
        q = "q{}".format(rid)
        lines = ["  const int {q} = rv{r} ? {pos} + ({off}) : {pos};".format(q=q, r=rid, pos=pos, off=off)]
        if lay.outer == "i" and dj:
            lines.append("  const int c{r} = rv{r} ? j + ({dj}) : j;".format(r=rid, dj=dj))
            rest = " + c{} * {}".format(rid, NK)
        lines.append("  const {ft}* __restrict__ p{r} = sf_cl_map({s} + ({q} - ({q} / {P}) * {P}) * {pl}{rest}, {q} / {P});"
                     .format(q=q, r=rid, ft=ft, s=slot, P=lay.P, pl=lay.plane, rest=rest))
        return "\n".join(lines)

    def _address(self, field, prow, kk):
        if field in self.layout.slot and self.layout.outer == "k":
            return "sf_cl_at<{}, {}, {}>({}, {})".format(
                ctype_of(self.program.fields[field].data_type), self.layout.P, self.layout.C, prow, kk)
        return super()._address(field, prow, kk)

    def _element(self, field, prow, kk):
        if field in self.layout.slot and self.layout.outer == "k":
            return "*" + self._address(field, prow, kk)
        return super()._element(field, prow, kk)


def generate(program, layout, specialize=None):
    """(kernel name, source, launch args) of the cluster kernel of ``program``."""
    fields = program.fields
    lay = layout
    T = lay.threads
    NI, NJ, NK = program.shape3
    gfields = lay.inputs + [o for o in program.outputs]
    gname = {f: "g{}".format(n) for n, f in enumerate(gfields)}
    scalars = []
    gens = []
    for op in program.ops:
        gen = ClusterOpGen(op, program, lay, specialize)
        gens.append(gen)
        scalars += [s for s in gen.scalars if s not in scalars]
    sname = {s: "sc{}".format(n) for n, s in enumerate(scalars)}
    params = ["const {}* __restrict__ {}".format(ctype_of(fields[f].data_type), gname[f]) for f in lay.inputs]
    params += ["{}* __restrict__ {}".format(ctype_of(fields[f].data_type), gname[f]) for f in program.outputs]
    params += ["const {} {}".format(ctype_of(fields[s].data_type), sname[s]) for s in scalars]

    body = ["  extern __shared__ __align__(16) unsigned char sf_smem[];",
            "  const int lo = (int)sf_cluster_rank() * {};".format(lay.P),
            "  const int n_own = min({}, lo + {}) - lo;".format(lay.n, lay.P)]
    sm = {f: "sm{}".format(n) for n, f in enumerate(lay.smem)}
    for f in lay.smem:
        ft = ctype_of(fields[f].data_type)
        body.append("  {}* const {} = reinterpret_cast<{}*>(sf_smem + {});".format(ft, sm[f], ft, lay.offset[f]))
    # full-dimensional inputs -> the owner's shared memory, 16-byte vectors where every range allows them
    for f in lay.loaded:
        ft, nb = ctype_of(fields[f].data_type), fields[f].data_type.bytes
        vl = max(1, 16 // nb)
        if (lay.P * lay.plane) % vl or (lay.n * lay.plane) % vl:
            vl = 1
        body.append("  for (int e = threadIdx.x * {vl}; e < n_own * {pl}; e += {step})\n"
                    "    *reinterpret_cast<SfVec<{ft}, {vl}>*>({s} + e) = "
                    "*reinterpret_cast<const SfVec<{ft}, {vl}>*>({g} + (i64)lo * {pl} + e);".format(
                        vl=vl, pl=lay.plane, step=T * vl, ft=ft, s=sm[f], g=gname[f]))
    for m, (op, gen) in enumerate(zip(program.ops, gens)):
        if m in lay.barriers:
            body.append("  sf_cluster_sync();")
        V = gen.V
        kv = NK // V
        body.append("  {{   // {}".format(op.name))
        for f in gen.in_fields:
            if f in gname and f not in lay.slot:
                body.append("  const {}* __restrict__ {} = {};".format(
                    ctype_of(fields[f].data_type), gen.canon[f], gname[f]))
        if op.name in gname:
            body.append("  {}* __restrict__ fout = {};".format(ctype_of(op.data_type), gname[op.name]))
        body.append("  for (int it = threadIdx.x; it < n_own * {} / {}; it += {}) {{".format(lay.plane, V, T))
        if lay.outer == "i":
            body.append("  const int k0 = (it % {}) * {}; const int j = (it / {}) % {}; const int i = lo + it / {};".format(
                kv, V, kv, NJ, kv * NJ))
        elif lay.outer == "j":
            body.append("  const int k0 = (it % {}) * {}; const int j = lo + it / {}; const int i = 0;".format(kv, V, kv))
        else:
            body.append("  const int k0 = lo + it * {}; const int j = 0; const int i = 0;".format(V))
        body.append("  (void)i; (void)j;")
        for s in gen.scalars:
            body.append("  const {} {} = sf_keep({});".format(ctype_of(fields[s].data_type), gen.scanon[s], sname[s]))
        cell, lines, results = gen.emit_cell()
        body += cell + lines + [gen.result_line(results)]
        ot = ctype_of(op.data_type)
        if op.name in lay.slot:
            body.append("  sf_stv<{}, {}>({} + it * {}, res);".format(ot, V, sm[op.name], V))
        if op.name in gname:
            body.append("  sf_stv<{}, {}>(fout + ({}), res);".format(ot, V, gen.out_index()))
        body.append("  }")
        body.append("  }")
    body.append("  sf_cluster_sync();          // no CTA leaves while a peer may still read its shared memory")
    text = "\n".join(body)
    digest = hashlib.sha1((text + ";".join(params) + repr((lay.C, T))).encode()).hexdigest()[:12]
    name = "sf_cluster_{}".format(digest)
    src = ('extern "C" __global__ void __cluster_dims__({}, 1, 1) __launch_bounds__({})\n{}({})\n{{\n{}\n}}\n'.format(
        lay.C, T, name, ", ".join(params), text))
    args = [("buf", f) for f in gfields] + [("scalar", fields[s].data_type, s) for s in scalars]
    return name, src, args


def lower_program_cluster(lowered, layout, specialize=None) -> LaunchSpec:
    """The whole program as one launch of one cluster (``layout.fits`` must hold)."""
    program = lowered.program
    name, src, args = generate(program, layout, specialize)
    block = (layout.threads, 1, 1)
    lowered.kernels[name] = KernelSpec(name, src, block, "cluster")
    C = layout.C
    launch = LaunchSpec(kernel=name, grid_fn=lambda b, e: (C, 1, 1), block=block, smem=layout.smem_bytes,
                        args=args, ops=[op.name for op in program.ops], reads=list(layout.inputs),
                        writes=list(program.outputs), cells_per_unit=program.cells, family="cluster",
                        info=layout.describe())
    lowered.launches.append(launch)
    return launch
